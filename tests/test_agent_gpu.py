"""End-to-end GPU parity: the B200 A2CAgent (CUDA kernels through the C ABI) vs
 (a) the committed golden fixtures produced by the REAL reference A2CAgent (tests/golden/agent_*.pt) and
 (b) the CPU oracle at a larger shape,
on identical env tapes, initial weights and sampling noise.  fp32 path (mixed_precision: False).

Tolerances: rollout tensors / normalised batch: rtol 1e-4; per-minibatch losses / KL: rtol 2e-3;
weights after 2 epochs (8-16 Adam steps): atol 2e-5 (Adam divides by sqrt(v): tiny-gradient elements
amplify 1e-7 differences); lr sequence and running-stat counts: exact.
"""
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as O

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')
DEV = 'cuda:0'
RUNS = tempfile.TemporaryDirectory(prefix='b200_test_runs_')      # the agents' train_dir: private to this process, removed at exit


class TapeEnvGPU:
    """GPU twin of oracle.ppo_oracle.TapeEnv / tests/golden/gen_golden.py::TapeVecEnv."""

    def __init__(self, obs_tape, done_tape, timeout_tape, A, autoreset='same_step', act_bounds=(-1.0, 1.0)):
        self.obs_tape, self.done_tape, self.timeout_tape = obs_tape.to(DEV), done_tape.to(DEV), timeout_tape.to(DEV)
        self.A, self.autoreset, self.i, self.act_bounds = A, autoreset, 0, act_bounds

    def reset(self):
        self.i = 0
        return self.obs_tape[0].clone()

    def step(self, actions):
        rew = -(actions * actions).sum(-1) * 0.1
        self.i += 1
        j = self.i % self.obs_tape.shape[0]
        return self.obs_tape[j].clone(), rew, self.done_tape[j].clone(), {'time_outs': self.timeout_tape[j].clone()}

    def get_env_info(self):
        from rl_games_b200.common import Box
        info = {'observation_space': Box(-np.inf, np.inf, (self.obs_tape.shape[-1],)), 'action_space': Box(self.act_bounds[0], self.act_bounds[1], (self.A,))}
        if self.autoreset != 'same_step':
            info['autoreset_mode'] = self.autoreset
        return info

    def get_env_state(self):
        return None

    def set_env_state(self, s):
        pass


def make_agent(cfg_over, N, H, D, A, units, mb, env, init_state, rnn_units=0, rnn_before_mlp=True, activation='elu', space_over=None, network_over=None):
    from rl_games_b200.runner import Runner
    network = {'name': 'actor_critic', 'separate': False,
               'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None', 'mu_init': {'name': 'default'},
                                        'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
               'mlp': {'units': list(units), 'activation': activation, 'initializer': {'name': 'default'}}}
    network['space']['continuous'].update(space_over or {})          # e.g. min_sigma (agent_minsigma.pt)
    network.update(network_over or {})                               # e.g. separate: True (agent_separate.pt)
    if rnn_units:
        network['rnn'] = {'name': 'lstm', 'units': rnn_units, 'layers': 1, 'before_mlp': rnn_before_mlp}
    config = {'name': 'gpu_parity', 'env_name': 'unused', 'reward_shaper': {'scale_value': 1.0}, 'device': DEV,
              'multi_gpu': False, 'mixed_precision': False, 'normalize_input': True, 'normalize_value': True,
              'value_bootstrap': True, 'normalize_advantage': True, 'gamma': 0.99, 'tau': 0.95, 'learning_rate': 3e-4,
              'lr_schedule': 'adaptive', 'kl_threshold': 0.008, 'grad_norm': 1.0, 'entropy_coef': 0.0, 'truncate_grads': True,
              'e_clip': 0.2, 'clip_value': True, 'use_smooth_clamp': True, 'bound_loss_type': 'regularisation',
              'bounds_loss_coef': 0.0, 'max_epochs': 100, 'num_actors': N, 'horizon_length': H, 'minibatch_size': mb,
              'mini_epochs': 4, 'critic_coef': 2, 'print_stats': False, 'train_dir': RUNS.name}
    config.update(cfg_over)
    config['env_info'] = env.get_env_info()
    config['vec_env'] = env
    params = {'seed': 7, 'algo': {'name': 'a2c_continuous'}, 'model': {'name': 'continuous_a2c_logstd'}, 'network': network,
              'config': config}
    r = Runner()
    r.load({'params': params})
    r.params['config']['vec_env'] = env
    agent = r.algo_factory.create(r.algo_name, base_name='parity', params=r.params)
    agent.model.load_state_dict({k: v.to(DEV) for k, v in init_state.items()}, strict=False)
    agent.init_tensors()
    agent._repack()
    agent.obs = agent.env_reset()
    return agent


def _check_epoch(agent, ref_state, ref_ds, ref_losses, ref_lr, units, tight=True, lstm=False):
    fl = O.swap_and_flatten01
    torch.testing.assert_close(fl(agent.advs_n).cpu(), ref_ds['advantages'], rtol=2e-4, atol=2e-5)
    torch.testing.assert_close(fl(agent.returns_n.unsqueeze(2)).cpu(), ref_ds['returns'], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(fl(agent.old_values_n.unsqueeze(2)).cpu(), ref_ds['old_values'], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(fl(agent.neglogpacs).cpu(), ref_ds['old_logp_actions'], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(fl(agent.actions).cpu(), ref_ds['actions'], rtol=1e-5, atol=1e-5)
    if ref_ds.get('rnn_masks') is not None:
        assert torch.equal(fl(agent.valid).cpu(), ref_ds['rnn_masks'])
    st = agent.last_stats
    for col, key in ((0, 'a'), (1, 'c'), (2, 'e'), (4, 'kl')):
        if ref_losses.get(key) is not None:
            torch.testing.assert_close(st[:, col], ref_losses[key], rtol=2e-3, atol=2e-6, msg=lambda m: key + ': ' + m)
    assert agent.last_lr == pytest.approx(ref_lr, rel=1e-12)
    sd = agent.model.state_dict()
    for k in O.param_names(len(units), lstm=lstm, separate=getattr(agent.model, 'separate', False)):
        torch.testing.assert_close(sd[k].cpu(), ref_state[k], rtol=1e-3, atol=2e-5, msg=lambda m: k + ': ' + m)
    for pre in ('running_mean_std.', 'value_mean_std.'):
        if pre + 'count' not in ref_state:          # that normaliser is switched off in this fixture: same key set as the reference
            assert pre + 'count' not in sd
            continue
        assert int(sd[pre + 'count']) == int(ref_state[pre + 'count'])
        torch.testing.assert_close(sd[pre + 'running_mean'].cpu(), ref_state[pre + 'running_mean'].reshape(-1), rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(sd[pre + 'running_var'].cpu(), ref_state[pre + 'running_var'].reshape(-1), rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize('name', ['agent_base.pt', 'agent_masked.pt', 'agent_hardclip.pt', 'agent_lstm.pt', 'agent_rmsadv.pt'])
@pytest.mark.parametrize('graph', [False, True])
def test_agent_matches_reference_golden(name, graph):
    _golden_run(name, graph)


@pytest.mark.parametrize('graph', [False, True])
def test_lstm_after_mlp_agent_matches_reference_golden(graph):
    """rnn before_mlp: False, the reference default (network_builder.py:253-272): same kernels as agent_lstm.pt, composed
    trunk -> LSTM window -> heads; the fixture comes from the reference itself (tests/golden/gen_golden.py lstm_after)"""
    _golden_run('agent_lstm_after.pt', graph, {})


@pytest.mark.parametrize('graph', [False, True])
def test_standard_schedule_agent_matches_reference_golden(graph):
    """schedule_type 'standard' (what the shipped mjlab configs use): the adaptive-KL scheduler steps once per mini-epoch on the mean
    KL, inside the optimiser kernel of the mini-epoch's last minibatch -- also when the update phase replays as a CUDA graph"""
    _golden_run('agent_sched_standard.pt', graph, {})


@pytest.mark.parametrize('name', ['agent_misc.pt', 'agent_rescale.pt', 'agent_minsigma.pt'])
@pytest.mark.parametrize('graph', [False, True])
def test_agent_matches_reference_golden_more_config_keys(name, graph):
    """agent_misc.pt: linear LR + entropy schedule (first minibatch of an epoch on the previous epoch's value), all normalisers off,
    full reward shaper, unclipped actions into a non-unit box; agent_rescale.pt: ppo: False, clip + rescale into that box, masked
    rows, bound loss; agent_minsigma.pt: the sigma floor of the 'exp' parametrisation (models.py:296-300; configs/mjlab/ppo_lift_cube_yam.yaml):
    the kernels read log(exp(raw) + min_sigma) and their log-std gradient is chained to the raw parameter, with an entropy bonus (whose
    gradient reaches only sigma), hard clip, bound loss, unclipped actions, masked rows.  Validated kernels, flag combinations no other
    GPU test sets."""
    _golden_run(name, graph)


@pytest.mark.parametrize('name', ['agent_lstm_masked.pt', 'agent_lstm_after_masked.pt'])
@pytest.mark.parametrize('graph', [False, True])
def test_lstm_on_next_step_autoreset_env_matches_reference_golden(name, graph):
    """envpool-style envs with an LSTM policy (a2c_common.py:1097-1106, :1180-1191): masked filler rows, the absorbed state re-zeroed in
    the rollout, the train-time reset also entering the first real row"""
    _golden_run(name, graph, {})


def _golden_run(name, graph, extra=None):
    g = torch.load(os.path.join(GOLDEN, name), weights_only=False)
    cfgk = g['config']
    over = {k: cfgk[k] for k in ('clip_value', 'use_smooth_clamp', 'bound_loss_type', 'bounds_loss_coef', 'entropy_coef',
                                 'truncate_grads', 'value_bootstrap', 'mini_epochs', 'lr_schedule', 'weight_decay', 'critic_coef', 'seq_length',
                                 'normalize_rms_advantage', 'adv_rms_momentum', 'schedule_type', 'learning_rate', 'kl_threshold',
                                 'max_epochs', 'schedule_entropy', 'normalize_input', 'normalize_value', 'normalize_advantage', 'clip_actions',
                                 'games_to_track', 'e_clip', 'tau', 'gamma', 'ppo')
            if k in cfgk}
    over.setdefault('lr_schedule', None)
    over['b200_cuda_graph'] = graph
    if g.get('reward_shaper'):
        over['reward_shaper'] = dict(g['reward_shaper'])
    over.update(extra or {})
    env = TapeEnvGPU(g['obs_tape'], g['done_tape'], g['timeout_tape'], g['A'], g['autoreset'], g.get('act_bounds', (-1.0, 1.0)))
    lstm = g.get('rnn_units', 0) > 0
    agent = make_agent(over, g['N'], g['H'], g['D'], g['A'], g['units'], g['mb'], env, g['init_state'], rnn_units=g.get('rnn_units', 0),
                       rnn_before_mlp=bool(g.get('rnn_before_mlp', True)), space_over=g.get('space_over'), network_over=g.get('network_over'))
    for ep, ref in enumerate(g['epochs_out']):
        agent.epoch_num += 1
        agent.train_epoch(noise=g['noise'][ep].to(DEV))
        assert torch.equal(agent.dones_buf.cpu(), ref['mb_dones'])
        torch.testing.assert_close(agent.rewards.cpu().unsqueeze(2), ref['mb_rewards'], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(agent.values.cpu().unsqueeze(2), ref['mb_values'], rtol=1e-4, atol=1e-5)
        nmb = agent.num_minibatches
        # reference returns per-minibatch a/c/entropy lists, per-mini-epoch mean KLs
        st = agent.last_stats
        torch.testing.assert_close(torch.stack([st[e * nmb:(e + 1) * nmb, 4].mean() for e in range(agent.mini_epochs_num)]),
                                   ref['kls'], rtol=2e-3, atol=2e-6)
        _check_epoch(agent, ref['state'], ref['dataset'], {'a': ref['a_losses'], 'c': ref['c_losses'], 'e': ref['entropies']},
                     ref['last_lr'], g['units'], lstm=lstm)
        torch.testing.assert_close(agent.game_rewards.mean, ref['game_rewards_mean'].reshape(-1), rtol=1e-4, atol=1e-5)
        assert agent.game_rewards.current_size == ref['game_rewards_size']
        torch.testing.assert_close(agent.game_lengths.mean, ref['game_lengths_mean'].reshape(-1), rtol=1e-5, atol=1e-5)
    return agent


@pytest.mark.parametrize('masked', [False, True])
def test_agent_matches_oracle_medium(masked):
    """N=256, H=16, D=60, A=8, MLP[64,32,16], mb=1024: exercises multi-block kernels and chunked minibatch rows."""
    N, H, D, A, units, mb, epochs = 256, 16, 60, 8, [64, 32, 16], 1024, 2
    obs_tape, done_tape, tout_tape = O.make_tapes(H * epochs + 1, N, D, seed=11)
    params = O.init_params(D, units, A, seed=3)
    g = torch.Generator().manual_seed(5)
    for k in params:
        if k.endswith('bias') or k.endswith('sigma'):
            params[k] = params[k] + torch.randn(params[k].shape, generator=g) * 0.05
    noise = torch.randn(epochs, H, N, A, generator=g)
    cfg = {'mask_autoreset_rows': masked, 'mini_epochs': 2}
    oag = O.OracleAgent(O.TapeEnv(obs_tape, done_tape, tout_tape), params, D, A, units, N, H, mb, cfg)
    oag.obs = oag.env_reset()
    env = TapeEnvGPU(obs_tape, done_tape, tout_tape, A, 'next_step' if masked else 'same_step')
    agent = make_agent({'mini_epochs': 2}, N, H, D, A, units, mb, env, params)
    for ep in range(epochs):
        out = oag.train_epoch(noise[ep])
        agent.epoch_num += 1
        agent.train_epoch(noise=noise[ep].to(DEV))
        ref_state = {k: v.detach() for k, v in oag.model.p.items()}
        for pre, m in (('running_mean_std.', oag.model.running_mean_std), ('value_mean_std.', oag.model.value_mean_std)):
            ref_state[pre + 'running_mean'], ref_state[pre + 'running_var'], ref_state[pre + 'count'] = \
                m.running_mean, m.running_var, m.count
        ds = {k: oag.dataset[k] for k in ('advantages', 'returns', 'old_values', 'old_logp_actions', 'actions', 'rnn_masks')}
        _check_epoch(agent, ref_state, ds, {'a': torch.stack(out['a_loss']), 'c': torch.stack(out['c_loss']),
                                            'e': torch.stack(out['entropy']), 'kl': torch.stack(out['kl'])}, oag.last_lr, units)


def test_checkpoint_roundtrip_and_reference_keys(tmp_path):
    N, H, D, A, units, mb = 64, 8, 6, 3, [16, 8], 128
    obs_tape, done_tape, tout_tape = O.make_tapes(H * 3 + 1, N, D, seed=2)
    env = TapeEnvGPU(obs_tape, done_tape, tout_tape, A)
    agent = make_agent({}, N, H, D, A, units, mb, env, O.init_params(D, units, A, seed=1))
    agent.epoch_num += 1
    agent.train_epoch()
    fn = str(tmp_path / 'ckpt')
    agent.save(fn)
    ck = torch.load(fn + '.pth', weights_only=False)
    # reference checkpoint layout: a2c_common.py:825-850 + state-dict keys (SURVEY 8b)
    assert set(['model', 'epoch', 'frame', 'optimizer', 'last_mean_rewards']).issubset(ck.keys())
    exp = set(O.param_names(len(units))) | {p + s for p in ('running_mean_std.', 'value_mean_std.')
                                             for s in ('running_mean', 'running_var', 'count')}
    assert set(ck['model'].keys()) == exp
    assert ck['model']['running_mean_std.count'].shape == () and ck['model']['running_mean_std.count'].dtype == torch.int64
    assert len(ck['optimizer']['state']) == 1 + 2 * len(units) + 4
    env2 = TapeEnvGPU(obs_tape, done_tape, tout_tape, A)
    agent2 = make_agent({}, N, H, D, A, units, mb, env2, O.init_params(D, units, A, seed=9))
    agent2.restore(fn + '.pth')
    assert torch.equal(agent2.model.flat, agent.model.flat)
    assert torch.equal(agent2.model.exp_avg, agent.model.exp_avg)
    # reference semantics (a2c_common.py:852-866): the optimizer comes back with its lr (held for the first step after the restore),
    # the agent's own last_lr is not part of a checkpoint
    assert agent2._resume_opt_lr == agent.last_lr and agent2.last_lr == 3e-4 and agent2.epoch_num == agent.epoch_num
    assert agent2.get_full_state_weights()['optimizer']['param_groups'][0]['lr'] == agent.last_lr
    torch.testing.assert_close(agent2.opt_state[1:4], agent.opt_state[1:4], rtol=1e-12, atol=0)      # step, beta1^step, beta2^step


def test_resume_from_a_reference_checkpoint_continues_like_the_reference():
    """tests/golden/gen_golden.py resume: a checkpoint of the REAL reference loaded into a fresh trainer, one more epoch -> where the
    reference's own fresh agent landed (weights, adaptive LR, Adam step count, normaliser statistics, epoch / frame)"""
    g = torch.load(os.path.join(GOLDEN, 'agent_resume.pt'), weights_only=False)
    ref, ck = g['resumed_epoch'], g['checkpoint']
    env = TapeEnvGPU(g['obs_tape'], g['done_tape'], g['timeout_tape'], g['A'])
    agent = make_agent({'weight_decay': g['config']['weight_decay'], 'lr_schedule': 'adaptive'}, g['N'], g['H'], g['D'], g['A'], g['units'], g['mb'],
                       env, g['init_state'])
    agent.set_full_state_weights({k: ({kk: vv.to(DEV) for kk, vv in v.items()} if k == 'model' else v) for k, v in ck.items()})
    agent.obs = agent.env_reset()
    agent.epoch_num += 1
    agent.train_epoch(noise=g['noise'][1].to(DEV))
    assert agent.epoch_num == ref['epoch_num'] and agent.frame == ref['frame']
    assert agent.last_lr == pytest.approx(ref['last_lr'], rel=1e-12)
    sd = agent.model.state_dict()
    for k in O.param_names(len(g['units'])):
        torch.testing.assert_close(sd[k].cpu(), ref['state'][k], rtol=1e-3, atol=2e-5, msg=lambda m: k + ': ' + m)
    out = agent.get_full_state_weights()
    assert float(out['optimizer']['state'][0]['step']) == ref['adam_step']


@pytest.mark.parametrize('mp', [False, True])
def test_masked_rows_contribute_zero_gradient(mp):
    """The reference's poison test (tests/test_ppo_masking.py:153-175), same call sequence: poison returns / values of the filler reset
    rows before prepare_dataset; one epoch of train_actor_critic from identical weights must give BIT-identical parameters (atol = 0) --
    masked value-normaliser moments, masked advantage normalisation, zero loss weight.  fp32 kernels and the bf16 tcgen05 kernels."""
    N, H, D, A, units, mb = (512, 8, 60, 8, [256, 128, 64], 2048) if mp else (64, 8, 6, 3, [16, 8], 128)
    obs_tape, done_tape, tout_tape = O.make_tapes(H + 1, N, D, seed=31)
    params = O.init_params(D, units, A, seed=5)
    g = torch.Generator().manual_seed(8)
    noise = torch.randn(H, N, A, generator=g).to(DEV)
    results = []
    for poison in (False, True):
        env = TapeEnvGPU(obs_tape, done_tape, tout_tape, A, autoreset='next_step')
        agent = make_agent({'mixed_precision': mp, 'mini_epochs': 2, 'b200_cuda_graph': False}, N, H, D, A, units, mb, env, params)
        # a first rollout so that the second one starts with pending reset rows at step 0 as well
        agent.play_steps(noise=noise)
        batch = agent.play_steps(noise=noise)
        garbage = batch['rnn_masks'] == 0.0
        assert 0 < int(garbage.sum()) < garbage.numel()
        if poison:
            batch['returns'] = batch['returns'].clone()
            batch['values'] = batch['values'].clone()
            batch['returns'][garbage] = 1e6
            batch['values'][garbage] = -1e6
        agent.set_train()
        agent.prepare_dataset(batch)
        for _ in range(agent.mini_epochs_num):
            for i in range(len(agent.dataset)):
                agent.train_actor_critic(agent.dataset[i])
        torch.cuda.synchronize()
        results.append({k: v.clone() for k, v in agent.model.state_dict().items()})
    clean, poisoned = results
    for k in clean:
        assert torch.equal(clean[k], poisoned[k]), f'parameter {k} differs: poisoned garbage rows leaked into the update'


def test_synthetic_env_training_runs_and_graph_replay_is_consistent():
    """c2-shaped (scaled down) synthetic env through the public Runner API; CUDA-graph replay vs eager updates
    from identical state must give identical weights (same kernels, same order => deterministic)."""
    from rl_games_b200.runner import Runner

    def build(graph):
        params = {'seed': 5, 'algo': {'name': 'a2c_continuous'}, 'model': {'name': 'continuous_a2c_logstd'},
                  'network': {'name': 'actor_critic', 'separate': False,
                              'space': {'continuous': {'mu_activation': 'None', 'sigma_activation': 'None',
                                                       'mu_init': {'name': 'default'},
                                                       'sigma_init': {'name': 'const_initializer', 'val': 0}, 'fixed_sigma': True}},
                              'mlp': {'units': [64, 32], 'activation': 'elu', 'initializer': {'name': 'default'}}},
                  'config': {'name': 'synt', 'env_name': 'b200_synthetic', 'reward_shaper': {'scale_value': 1.0}, 'device': DEV,
                             'normalize_input': True, 'normalize_value': True, 'normalize_advantage': True, 'gamma': 0.99,
                             'tau': 0.95, 'learning_rate': 3e-4, 'lr_schedule': 'adaptive', 'kl_threshold': 0.008,
                             'grad_norm': 1.0, 'entropy_coef': 0.0, 'truncate_grads': True, 'e_clip': 0.2, 'clip_value': True,
                             'use_smooth_clamp': True, 'bound_loss_type': 'regularisation', 'bounds_loss_coef': 0.0,
                             'num_actors': 1024, 'horizon_length': 16, 'minibatch_size': 4096, 'mini_epochs': 2,
                             'critic_coef': 2, 'print_stats': False, 'train_dir': RUNS.name,
                             'mixed_precision': False, 'b200_cuda_graph': graph,
                             'env_config': {'obs_dim': 60, 'act_dim': 8, 'device': DEV}}}
        r = Runner()
        r.load({'params': params})
        a = r.algo_factory.create(r.algo_name, base_name='synt', params=r.params)
        a.init_tensors()
        a.obs = a.env_reset()
        return a
    a, b = build(True), build(False)
    b.model.load_state_dict(a.model.state_dict())
    for _ in range(4):
        a.epoch_num += 1; b.epoch_num += 1
        a.train_epoch(); b.train_epoch()
    assert (a._graph_epoch is not None or a._graph_update is not None) and b._graph_update is None and b._graph_epoch is None
    assert torch.equal(a.model.flat, b.model.flat)
    assert a.last_lr == b.last_lr
    assert torch.isfinite(a.model.flat).all()
    assert a.game_rewards.current_size > 0


def test_bf16_tcgen05_agent_tracks_fp32_agent():
    """mixed_precision: True (bf16 tcgen05 kernels) vs mixed_precision: False (fp32 kernels) on the c2 architecture
    (obs 60, MLP [256,128,64], 8 actions), same tapes / weights / noise.  bf16 tolerance class (8-bit mantissa operands,
    fp32 accumulate): rollout outputs atol 5e-2, per-minibatch losses rtol 0.1 (+ small atol), parameter update
    direction cosine > 0.8 after one epoch of Adam steps."""
    _bf16_vs_fp32_agents(60, {})


@pytest.mark.parametrize('D', [256, 105])
def test_bf16_tcgen05_wide_agent_tracks_fp32_agent(D):
    """the same comparison on BASELINE configs[4]'s observation width (256) and a ragged one: layer 1 in its own kernels"""
    _bf16_vs_fp32_agents(D, {})


@pytest.mark.parametrize('extra', [{'ppo': False}, {'normalize_input': False, 'normalize_value': False, 'normalize_advantage': False},
                                   {'clip_actions': False}, {'clip_value': False, 'use_smooth_clamp': False},
                                   {'bounds_loss_coef': 0.001, 'bound_loss_type': 'bound'}, {'bounds_loss_coef': None},
                                   {'truncate_grads': False, 'weight_decay': 0.01, 'entropy_coef': 0.01}],
                         ids=lambda e: ','.join(f'{k}={v}' for k, v in e.items()))
def test_bf16_tcgen05_agent_tracks_fp32_agent_flag_matrix(extra):
    """every loss / shaping / optimiser flag the fused tcgen05 kernels branch on, against the fp32 kernels (which the reference golden
    runs pin): same tolerance class as the default comparison"""
    _bf16_vs_fp32_agents(60, dict(extra))


@pytest.mark.parametrize('D,units,activation', [(17, [128, 64, 32], 'relu'), (60, [128, 64, 32], 'tanh'), (111, [200, 100, 50], 'elu'), (60, [256, 128, 64], 'relu')])
def test_bf16_tcgen05_agent_other_geometries_and_activations_track_fp32_agent(D, units, activation):
    """three-layer MLPs narrower than the compiled tiles (zero-padded; [128, 64, 32] is configs/mujoco/walker2d.yaml) and relu / tanh
    networks on the tcgen05 kernels vs the fp32 kernels: the same tolerance class as the native geometry"""
    _bf16_vs_fp32_agents(D, {}, units=units, activation=activation)


def _bf16_vs_fp32_agents(D, extra, units=(256, 128, 64), activation='elu'):
    N, H, A, mb = 512, 8, 8, 2048
    units = list(units)
    obs_tape, done_tape, tout_tape = O.make_tapes(H + 1, N, D, seed=21)
    params = O.init_params(D, units, A, seed=4)
    g = torch.Generator().manual_seed(6)
    noise = torch.randn(H, N, A, generator=g).to(DEV)
    agents = []
    for mp in (False, True):
        env = TapeEnvGPU(obs_tape, done_tape, tout_tape, A)
        a = make_agent({'mixed_precision': mp, 'mini_epochs': 2, 'b200_cuda_graph': False, **extra}, N, H, D, A, units, mb, env, params, activation=activation)
        assert a.use_tc == mp and getattr(a, 'tc_wide', False) == (mp and D > 64)
        a.epoch_num += 1
        a.train_epoch(noise=noise)
        agents.append(a)
    f, t = agents
    torch.testing.assert_close(t.values, f.values, rtol=0, atol=6e-2)
    torch.testing.assert_close(t.mus, f.mus, rtol=0, atol=6e-2)   # after the update: last mini-epoch's mu write-back
    torch.testing.assert_close(t.advs_n, f.advs_n, rtol=0, atol=0.15)
    sf, st = f.last_stats, t.last_stats
    torch.testing.assert_close(st[:, 0], sf[:, 0], rtol=0.1, atol=2e-2)     # a_loss
    torch.testing.assert_close(st[:, 1], sf[:, 1], rtol=0.1, atol=2e-2)     # c_loss
    torch.testing.assert_close(st[:, 2], sf[:, 2], rtol=1e-3, atol=1e-3)    # entropy (depends on sigma only)
    torch.testing.assert_close(st[:, 4], sf[:, 4], rtol=0.35, atol=3e-4)    # kl
    init = torch.cat([params[k].reshape(-1) for k in O.param_names(3)])
    # flat order differs from param_names order only by the head packing; compare per tensor through state_dict
    sdf, sdt = f.model.state_dict(), t.model.state_dict()
    for k in O.param_names(3):
        if k.endswith('weight'):
            du_f = (sdf[k].cpu() - params[k]).flatten(); du_t = (sdt[k].cpu() - params[k]).flatten()
            cos = float(du_f @ du_t / (du_f.norm() * du_t.norm() + 1e-20))
            assert cos > 0.8, (k, cos)
    assert 0.4 < t.last_lr / f.last_lr < 2.5
    if t.normalize_input:
        assert int(t.model.running_mean_std.count) == int(f.model.running_mean_std.count)


@pytest.mark.parametrize('opt', [{'b200_pdl': True}, {'b200_pipelined_wgrad': True}, {'b200_pdl': True, 'b200_cuda_graph': True}])
def test_tc_agent_launch_options_do_not_change_results(opt):
    """programmatic dependent launch (b200_pdl) only changes WHEN the chain kernels may start, never what they compute: weights
    after two epochs are bit-identical to the plain stream-ordered run (eager and whole-epoch graph).  The pipelined
    weight-gradient kernel (b200_pipelined_wgrad) sums rows in 64-row halves: fp32 accumulation-order agreement."""
    from rl_games_b200 import ops
    N, H, D, A, units, mb = 1024, 8, 60, 8, [256, 128, 64], 4096
    obs_tape, done_tape, tout_tape = O.make_tapes(2 * H + 1, N, D, seed=23)
    params = O.init_params(D, units, A, seed=5)
    g = torch.Generator().manual_seed(7)
    noise = [torch.randn(H, N, A, generator=g).to(DEV) for _ in range(2)]
    out = []
    try:
        for over in ({}, opt):
            env = TapeEnvGPU(obs_tape, done_tape, tout_tape, A)
            cfg = {'mixed_precision': True, 'mini_epochs': 2, 'b200_cuda_graph': False}
            cfg.update(over)
            a = make_agent(cfg, N, H, D, A, units, mb, env, params)
            assert a.use_tc
            for e in range(2):
                a.epoch_num += 1
                a.train_epoch(noise=noise[e])
            torch.cuda.synchronize()
            out.append((a.model.flat.clone(), a.last_stats.clone(), a.last_lr))
    finally:
        ops.set_pdl(False)
    (f0, s0, lr0), (f1, s1, lr1) = out
    assert torch.isfinite(f1).all()
    if 'b200_pipelined_wgrad' in opt:
        torch.testing.assert_close(f1, f0, rtol=0, atol=2e-4)        # Adam steps of 3e-4: a sign flip of a ~0 gradient moves a weight by <= lr
        torch.testing.assert_close(s1[:, :5], s0[:, :5], rtol=2e-2, atol=1e-3)
    else:
        assert torch.equal(f1, f0) and torch.equal(s1, s0) and lr1 == lr0


@pytest.mark.parametrize('name,N,H,D,A,mb,masked,mp', [
    ('c3_ant_envpool_shape', 4096, 64, 27, 8, 32768, True, False),     # BASELINE configs[2]: next_step autoreset => masked path
    ('c5_per_gpu_shape', 16384, 32, 256, 8, 32768, False, False),      # BASELINE configs[4] per-GPU shard (obs 256): fp32 path
    ('c2_shape_bf16', 16384, 16, 60, 8, 32768, False, True),           # BASELINE configs[1] on the tcgen05 path
])
def test_full_size_configs_one_epoch_vs_oracle(name, N, H, D, A, mb, masked, mp):
    """BASELINE.json full-size shapes: one complete epoch (rollout -> GAE -> 1 mini-epoch of updates) against the CPU oracle
    on identical tapes / weights / noise.  fp32 path: rollout + normalised batch rtol 1e-4, losses rtol 5e-3, weights atol 5e-5;
    bf16 path: bf16 tolerance class."""
    units = [256, 128, 64]
    g = torch.Generator().manual_seed(17)
    T = H + 1
    obs_tape = torch.randn(T, N, D, generator=g) * 1.5 + 0.3
    done_tape = (torch.rand(T, N, generator=g) < 0.03).to(torch.uint8)
    tout_tape = (torch.rand(T, N, generator=g) < 0.3) & done_tape.bool()
    params = O.init_params(D, units, A, seed=6)
    noise = torch.randn(H, N, A, generator=g)
    oag = O.OracleAgent(O.TapeEnv(obs_tape, done_tape, tout_tape), params, D, A, units, N, H, mb,
                        {'mask_autoreset_rows': masked, 'mini_epochs': 1}, matmul_dtype=torch.bfloat16 if mp else None)
    oag.obs = oag.env_reset()
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    out = oag.train_epoch(noise)
    env = TapeEnvGPU(obs_tape, done_tape, tout_tape, A, 'next_step' if masked else 'same_step')
    agent = make_agent({'mini_epochs': 1, 'mixed_precision': mp}, N, H, D, A, units, mb, env, params)
    agent.epoch_num += 1
    agent.train_epoch(noise=noise.to(DEV))
    fl = O.swap_and_flatten01
    st = agent.last_stats
    if not mp:
        assert torch.equal(agent.dones_buf.cpu(), oag.buf['dones'])
        torch.testing.assert_close(agent.values.cpu(), oag.buf['values'].squeeze(2), rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(fl(agent.advs_n).cpu(), oag.dataset['advantages'], rtol=1e-3, atol=1e-4)
        torch.testing.assert_close(st[:, 0], torch.stack(out['a_loss']), rtol=5e-3, atol=1e-5)
        torch.testing.assert_close(st[:, 1], torch.stack(out['c_loss']), rtol=5e-3, atol=1e-5)
        torch.testing.assert_close(st[:, 4], torch.stack(out['kl']), rtol=1e-2, atol=1e-6)
        assert agent.last_lr == pytest.approx(oag.last_lr, rel=1e-12)
        sd = agent.model.state_dict()
        for k in O.param_names(3):
            torch.testing.assert_close(sd[k].cpu(), oag.model.p[k].detach(), rtol=1e-3, atol=5e-5, msg=lambda m: k + ': ' + m)
        assert int(sd['running_mean_std.count']) == int(oag.model.running_mean_std.count)
        torch.testing.assert_close(sd['running_mean_std.running_mean'].cpu(), oag.model.running_mean_std.running_mean, rtol=1e-5, atol=1e-6)
    else:
        torch.testing.assert_close(agent.values.cpu(), oag.buf['values'].squeeze(2), rtol=0, atol=8e-2)
        torch.testing.assert_close(st[:, 0], torch.stack(out['a_loss']), rtol=0.15, atol=3e-3)
        torch.testing.assert_close(st[:, 1], torch.stack(out['c_loss']), rtol=0.1, atol=2e-2)
        torch.testing.assert_close(st[:, 4], torch.stack(out['kl']), rtol=0.3, atol=2e-4)
        assert int(agent.model.running_mean_std.count) == int(oag.model.running_mean_std.count)


def test_lstm_agent_matches_oracle_medium():
    """LSTM-before-MLP policy (BASELINE configs[3] structure, scaled down): N=128 envs, H=16, seq_length=4, obs 44, 5 actions, LSTM 32,
    MLP [64,32]; two epochs with episode ends inside the BPTT windows; fp32 path vs the CPU oracle (pinned to the reference by
    tests/golden/agent_lstm.pt)."""
    N, H, D, A, units, mb, hid, epochs = 128, 16, 44, 5, [64, 32], 512, 32, 2
    obs_tape, done_tape, tout_tape = O.make_tapes(H * epochs + 1, N, D, seed=31, p_done=0.08)
    params = O.init_params(D, units, A, seed=3, rnn_units=hid)
    g = torch.Generator().manual_seed(15)
    noise = torch.randn(epochs, H, N, A, generator=g)
    cfg = {'mini_epochs': 2, 'rnn_units': hid, 'seq_length': 4}
    oag = O.OracleAgent(O.TapeEnv(obs_tape, done_tape, tout_tape), params, D, A, units, N, H, mb, cfg)
    oag.obs = oag.env_reset()
    env = TapeEnvGPU(obs_tape, done_tape, tout_tape, A)
    agent = make_agent({'mini_epochs': 2, 'seq_length': 4}, N, H, D, A, units, mb, env, params, rnn_units=hid)
    assert agent.is_rnn and not agent.use_tc
    for ep in range(epochs):
        out = oag.train_epoch(noise[ep])
        agent.epoch_num += 1
        agent.train_epoch(noise=noise[ep].to(DEV))
        ref_state = {k: v.detach() for k, v in oag.model.p.items()}
        for pre, m in (('running_mean_std.', oag.model.running_mean_std), ('value_mean_std.', oag.model.value_mean_std)):
            ref_state[pre + 'running_mean'], ref_state[pre + 'running_var'], ref_state[pre + 'count'] = \
                m.running_mean, m.running_var, m.count
        ds = {k: oag.dataset[k] for k in ('advantages', 'returns', 'old_values', 'old_logp_actions', 'actions', 'rnn_masks')}
        _check_epoch(agent, ref_state, ds, {'a': torch.stack(out['a_loss']), 'c': torch.stack(out['c_loss']),
                                            'e': torch.stack(out['entropy']), 'kl': torch.stack(out['kl'])}, oag.last_lr, units, lstm=True)
        # rollout-side state snapshots (mb_rnn_states, a2c_common.py:1081-1083) and the carried states
        torch.testing.assert_close(agent.rnn_h0.cpu(), oag.mb_rnn_states[0].squeeze(1), rtol=1e-4, atol=1e-5)
        torch.testing.assert_close(agent.rnn_c0.cpu(), oag.mb_rnn_states[1].squeeze(1), rtol=1e-4, atol=1e-5)
        torch.testing.assert_close(agent.rnn_h.cpu(), oag.rnn_states[0][0], rtol=1e-4, atol=1e-5)


def test_lstm_c4_geometry_full_width_vs_oracle():
    """BASELINE configs[3] geometry at full width: 8192 envs, obs 348, 17 actions (Humanoid-v5), LSTM 256 before the MLP [512, 256, 128]
    (configs/mujoco/humanoid_envpool.yaml:23), seq_length 4 -- horizon 8 (two BPTT windows per env; the horizon only repeats windows), one
    mini-epoch of 4 minibatches, fp32 kernels vs the CPU oracle on identical tapes / weights / noise: rollout values and states rtol 1e-4,
    losses rtol 5e-3, weights atol 5e-5."""
    N, H, D, A, units, mb, hid = 8192, 8, 348, 17, [512, 256, 128], 16384, 256
    g = torch.Generator().manual_seed(41)
    T = H + 1
    obs_tape = torch.randn(T, N, D, generator=g) * 1.5 + 0.3
    done_tape = (torch.rand(T, N, generator=g) < 0.05).to(torch.uint8)
    tout_tape = (torch.rand(T, N, generator=g) < 0.3) & done_tape.bool()
    params = O.init_params(D, units, A, seed=9, rnn_units=hid)
    noise = torch.randn(H, N, A, generator=g)
    cfg = {'mini_epochs': 1, 'rnn_units': hid, 'seq_length': 4}
    oag = O.OracleAgent(O.TapeEnv(obs_tape, done_tape, tout_tape), params, D, A, units, N, H, mb, cfg)
    oag.obs = oag.env_reset()
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    out = oag.train_epoch(noise)
    env = TapeEnvGPU(obs_tape, done_tape, tout_tape, A)
    agent = make_agent({'mini_epochs': 1, 'seq_length': 4}, N, H, D, A, units, mb, env, params, rnn_units=hid)
    assert agent.is_rnn and not agent.use_tc and agent.model.rnn_units == hid
    agent.epoch_num += 1
    agent.train_epoch(noise=noise.to(DEV))
    st = agent.last_stats
    torch.testing.assert_close(agent.values.cpu(), oag.buf['values'].squeeze(2), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(agent.rnn_h.cpu(), oag.rnn_states[0][0], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(st[:, 0], torch.stack(out['a_loss']), rtol=5e-3, atol=1e-5)
    torch.testing.assert_close(st[:, 1], torch.stack(out['c_loss']), rtol=5e-3, atol=1e-5)
    torch.testing.assert_close(st[:, 4], torch.stack(out['kl']), rtol=1e-2, atol=1e-6)
    assert agent.last_lr == pytest.approx(oag.last_lr, rel=1e-12)
    sd = agent.model.state_dict()
    for k in O.param_names(3, lstm=True):
        torch.testing.assert_close(sd[k].cpu(), oag.model.p[k].detach(), rtol=1e-3, atol=5e-5, msg=lambda m: k + ': ' + m)


def test_rollout_precision_option_reproduces_the_fp32_rollout_exactly():
    """b200_rollout_fp32 (the reference's precision split: rollout outside autocast, a2c_common.py:581-600; update in bf16,
    a2c_continuous.py:173): with it the tcgen05 agent's rollout arena is BIT-identical to the fp32 agent's on the same weights / noise;
    without it (default: bf16 rollout, self-consistent with the bf16 update) the arena differs by the bf16 tolerance class, measured
    here: |dvalue| <= 6e-2, |dmu| <= 6e-2, and the first-minibatch importance ratio is exactly 1 only in the default mode."""
    N, H, D, A, units, mb = 512, 8, 60, 8, [256, 128, 64], 2048
    obs_tape, done_tape, tout_tape = O.make_tapes(H + 1, N, D, seed=33)
    params = O.init_params(D, units, A, seed=8)
    g = torch.Generator().manual_seed(9)
    noise = torch.randn(H, N, A, generator=g).to(DEV)
    ag = {}
    for name, cfg in (('fp32', {'mixed_precision': False}), ('tc', {'mixed_precision': True}),
                      ('tc_rollout_fp32', {'mixed_precision': True, 'b200_rollout_fp32': True})):
        # normalize_input off: the obs normaliser moves between the rollout and the first minibatch (model.train()), which would hide the precision effect
        a = make_agent({'mini_epochs': 1, 'b200_cuda_graph': False, 'normalize_input': False, **cfg}, N, H, D, A, units, mb,
                       TapeEnvGPU(obs_tape, done_tape, tout_tape, A), params)
        a._rollout(noise)
        a._gae_and_prepare()
        torch.cuda.synchronize()
        ag[name] = a
    f, t, tf = ag['fp32'], ag['tc'], ag['tc_rollout_fp32']
    assert tf.use_tc and tf.rollout_fp32 and not t.rollout_fp32
    for k in ('values', 'mus', 'neglogpacs', 'actions', 'rewards', 'advs_n', 'returns_n'):
        assert torch.equal(getattr(tf, k), getattr(f, k)), k
    torch.testing.assert_close(t.values, f.values, rtol=0, atol=6e-2)
    torch.testing.assert_close(t.mus, f.mus, rtol=0, atol=6e-2)
    # first minibatch: ratio = exp(old_neglogp - neglogp) == 1 <=> a_loss == -mean(adv) ... measured through the KL statistic (0 iff mu, sigma match)
    for a in (t, tf):
        a._minibatch_update(0, 0)
    torch.cuda.synchronize()
    kl_default, kl_split = float(t.stats[0, 4]), float(tf.stats[0, 4])
    # policy_kl of two IDENTICAL Gaussians is not 0 but A * (log(1 + 1e-5) + 1 / (2 (1 + 1e-5)) - 1/2) (the 1e-5 terms of torch_ext.py:27-36), sigma = 1 here
    import math
    kl_same = A * (math.log1p(1e-5) + 0.5 / (1.0 + 1e-5) - 0.5)
    assert abs(kl_default - kl_same) < 2e-6, (kl_default, kl_same)      # same arithmetic in rollout and update: the policy has not moved yet
    assert kl_default < kl_split < 5e-3, (kl_default, kl_split)          # fp32 behaviour policy vs bf16 re-evaluation: bf16 noise shows up as a spurious KL
    print('rollout precision: first-minibatch KL default (bf16 rollout) %.3e, reference split (fp32 rollout) %.3e' % (kl_default, kl_split))


@pytest.mark.parametrize('case', ['lstm_before_mlp', 'lstm_after_mlp', 'mlp_512_256_128', 'mlp_128_64_32_min_sigma'])
def test_layerwise_tensor_core_path_tracks_fp32_agent(case):
    """mixed_precision: True on an LSTM policy / an MLP wider than the fused tiles: every GEMM on the tensor cores (gemm_tc.cu, bf16
    operands, fp32 accumulate), the same host composition as the fp32 path.  Against the fp32 kernels on the same tapes / weights /
    noise: bf16 tolerance class (rollout outputs atol 6e-2, per-minibatch losses rtol 0.1, update direction cosine > 0.8).
    mlp_128_64_32_min_sigma: a geometry the FUSED kernels have, with a sigma floor (min_sigma; the fused kernels read the raw parameter from
    the packed arena, so the floored policy is routed layer by layer) -- the floor, its gradient chain and an entropy bonus on both paths."""
    N, H, D, A, mb = 256, 8, 44, 5, 1024
    units, rnn, before = ([64, 32], 32, True) if case == 'lstm_before_mlp' else (([64, 32], 32, False) if case == 'lstm_after_mlp' else ([512, 256, 128], 0, True))
    space_over, extra = None, {}
    if case == 'mlp_128_64_32_min_sigma':
        units, space_over, extra = [128, 64, 32], {'min_sigma': 0.2}, {'entropy_coef': 0.01}
    obs_tape, done_tape, tout_tape = O.make_tapes(H + 1, N, D, seed=51, p_done=0.08)
    params = O.init_params(D, units, A, seed=6, rnn_units=rnn, rnn_before_mlp=before)
    g = torch.Generator().manual_seed(16)
    noise = torch.randn(H, N, A, generator=g).to(DEV)
    agents = []
    for mp in (False, True):
        a = make_agent(dict({'mixed_precision': mp, 'mini_epochs': 2, 'b200_cuda_graph': False, 'seq_length': 4}, **extra), N, H, D, A, units, mb,
                       TapeEnvGPU(obs_tape, done_tape, tout_tape, A), params, rnn_units=rnn, rnn_before_mlp=before, space_over=space_over)
        assert a.gemm_tc == mp and not a.use_tc and a.model.min_sigma == (space_over or {}).get('min_sigma', 0.0)
        a.epoch_num += 1
        a.train_epoch(noise=noise)
        agents.append(a)
    f, t = agents
    torch.testing.assert_close(t.values, f.values, rtol=0, atol=6e-2)
    torch.testing.assert_close(t.mus, f.mus, rtol=0, atol=6e-2)
    sf, st = f.last_stats, t.last_stats
    torch.testing.assert_close(st[:, 0], sf[:, 0], rtol=0.1, atol=2e-2)
    torch.testing.assert_close(st[:, 1], sf[:, 1], rtol=0.1, atol=2e-2)
    torch.testing.assert_close(st[:, 4], sf[:, 4], rtol=0.35, atol=3e-4)
    sdf, sdt = f.model.state_dict(), t.model.state_dict()
    for k in O.param_names(len(units), lstm=bool(rnn)):
        if k.endswith('weight') or 'weight_' in k:
            du_f = (sdf[k].cpu() - params[k]).flatten(); du_t = (sdt[k].cpu() - params[k]).flatten()
            cos = float(du_f @ du_t / (du_f.norm() * du_t.norm() + 1e-20))
            assert cos > 0.8, (k, cos)
    if space_over:          # the floored sigma: the stored sigmas (rewritten by the last mini-epoch, datasets.py:33-43) are exp(raw) + min_sigma on
        # both paths -- equal up to what the two paths' slightly different updates did to raw (measured: 2e-6) -- and raw moved the same way
        torch.testing.assert_close(t.sigmas, f.sigmas, rtol=0, atol=1e-3)
        assert float(f.sigmas.min()) > space_over['min_sigma']
        ds_f, ds_t = sdf['a2c_network.sigma'].cpu() - params['a2c_network.sigma'], sdt['a2c_network.sigma'].cpu() - params['a2c_network.sigma']
        assert float(ds_f @ ds_t / (ds_f.norm() * ds_t.norm() + 1e-20)) > 0.8
